"""CUDA backend: drives the native sm_100a core for tensors that live on the GPU.

This is the layer the reference implements in mpi_xla_bridge_cuda.cpp (882 lines of
host C++ that synchronise the stream and hand pointers to MPI).  Here a communicator
owns peer-mapped HBM:

* a *control segment* (barrier flags, p2p rings, LL buffers, halo buffers) and
* a growable *staging segment* (+ its NVLS multicast alias),

both created with the CUDA VMM API inside ``libb2mpi.so``; the POSIX file descriptors
that name the physical allocations are exchanged between the local ranks over unix
domain sockets (``SCM_RIGHTS``), everything else over the gloo control plane.  Every
op is a kernel launch on the caller's current stream: nothing here synchronises the
host, so ops can be recorded into CUDA graphs (``mpi4jax_b200.jit``).
"""

from __future__ import annotations

import ctypes
import functools
import os
import socket
import sys
import tempfile
import threading
import uuid
import weakref
from typing import Optional

import torch
import torch.distributed as dist

from .. import native
from ..comm import ANY_SOURCE, ANY_TAG, Comm, MPIError, Status
from ..decorators import env_flag, env_float, env_int, setup_cuda_mpi
from ..native import codes

_MIN_STAGE = 64 << 20
_POISON = env_flag("MPI4JAX_B200_POISON", False)


class _RawDeviceBytes:
    """``__cuda_array_interface__`` view of raw device memory (for the poison debug mode)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False),
                                         "version": 2}


def _lib():
    if not native.HAS_CUDA_EXT:
        raise ImportError(
            "mpi4jax_b200: CUDA tensors need the native library, which failed to load "
            f"({native.CUDA_EXT_ERROR}); build it with `python -m mpi4jax_b200._src.native.build`."
        )
    return native.lib


def abort_or_raise(message: str, code: int = 1):
    """The reference's fail-fast path (mpi_ops_common.h:60-78): print
    ``r<rank> | MPI_<op> returned error code ... - aborting`` and kill the job."""
    sys.stderr.write(message + "\n")
    sys.stderr.flush()
    if env_flag("MPI4JAX_B200_ABORT_ON_ERROR", True):
        os._exit(code if 0 < code < 256 else 1)
    raise MPIError(message)


# ---------------------------------------------------------------------------
# control-plane helpers
# ---------------------------------------------------------------------------
def _all_gather_obj(comm: Comm, obj):
    out = [None] * comm.size
    if comm.size == 1:
        return [obj]
    dist.all_gather_object(out, obj, group=comm._group)
    return comm._in_rank_order(out)


def _exchange_fds(comm: Comm, fd: Optional[int]) -> dict:
    """Every rank that passes an fd sends a duplicate of it to all other ranks.
    Returns {source_rank: received_fd}."""
    if comm.size == 1:
        return {}
    token = uuid.uuid4().hex[:12]
    path = os.path.join(tempfile.gettempdir(), f"b2mpi-{os.getpid()}-{token}.sock")
    listener = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
    listener.bind(path)
    listener.listen(comm.size)
    info = _all_gather_obj(comm, (path, fd is not None))
    senders = [r for r, (_, has) in enumerate(info) if has and r != comm.rank]
    received: dict = {}
    errors: list = []

    def accept_all():
        try:
            for _ in senders:
                conn, _addr = listener.accept()
                with conn:
                    msg, fds, _flags, _a = socket.recv_fds(conn, 64, 1)
                    received[int(msg.decode())] = fds[0]
        except Exception as exc:  # pragma: no cover
            errors.append(exc)

    th = threading.Thread(target=accept_all, daemon=True)
    th.start()
    if fd is not None:
        for r, (peer_path, _) in enumerate(info):
            if r == comm.rank:
                continue
            with socket.socket(socket.AF_UNIX, socket.SOCK_STREAM) as s:
                s.connect(peer_path)
                socket.send_fds(s, [str(comm.rank).encode()], [fd])
    th.join(timeout=120)
    listener.close()
    try:
        os.unlink(path)
    except OSError:
        pass
    if errors or th.is_alive():
        raise MPIError(f"file-descriptor exchange failed: {errors}")
    dist.barrier(group=comm._group)
    return received


class _Segment:
    """A symmetric segment (+ optional multicast alias) shared by all ranks of a comm."""

    def __init__(self, comm: Comm, device: int, nbytes: int, mode: str, want_mc: bool):
        lib = _lib()
        self.comm = comm
        self.seg = None
        self.mc = None
        mode_code = 0 if mode == "vmm" else 1
        seg = lib.b2_seg_create(device, comm.rank, comm.size, nbytes, mode_code)
        oks = _all_gather_obj(comm, bool(seg))
        if not all(oks):
            err = native.last_error()
            if seg:
                lib.b2_seg_destroy(seg)
            raise MPIError(f"symmetric segment allocation failed on ranks "
                           f"{[r for r, ok in enumerate(oks) if not ok]}: {err}")
        self.seg = seg
        self.bytes = int(lib.b2_seg_bytes(seg))
        if comm.size > 1:
            if mode == "vmm":
                fd = lib.b2_seg_export_fd(seg)
                if fd < 0:
                    raise MPIError(f"exporting the segment failed: {native.last_error()}")
                for peer, pfd in _exchange_fds(comm, fd).items():
                    rc = lib.b2_seg_import_fd(seg, peer, pfd)
                    os.close(pfd)
                    if rc != 0:
                        raise MPIError(f"mapping rank {peer}'s segment failed: {native.last_error()}")
            else:
                buf = ctypes.create_string_buffer(64)
                if lib.b2_seg_ipc_handle(seg, buf) != 0:
                    raise MPIError(f"cudaIpcGetMemHandle failed: {native.last_error()}")
                handles = _all_gather_obj(comm, bytes(buf.raw))
                for peer, h in enumerate(handles):
                    if peer == comm.rank:
                        continue
                    hb = ctypes.create_string_buffer(h, 64)
                    if lib.b2_seg_import_ipc(seg, peer, hb) != 0:
                        raise MPIError(f"cudaIpcOpenMemHandle failed: {native.last_error()}")
            dist.barrier(group=comm._group)
        if want_mc and mode == "vmm" and comm.size > 1:
            self._setup_multicast(device)

    def _setup_multicast(self, device: int) -> None:
        lib = _lib()
        comm = self.comm
        mc = None
        fd = None
        if comm.rank == 0:
            mc = lib.b2_mc_create(device, comm.size, self.bytes)
            if mc:
                fd = lib.b2_mc_export_fd(mc)
                if fd < 0:
                    lib.b2_mc_destroy(mc)
                    mc, fd = None, None
        ok0 = _all_gather_obj(comm, bool(mc) if comm.rank == 0 else True)[0]
        if not ok0:
            return                      # multicast unavailable: plain P2P paths only
        got = _exchange_fds(comm, fd)
        if comm.rank != 0:
            mc = lib.b2_mc_import(device, got[0], self.bytes)
            os.close(got[0])
        ok = bool(mc) and lib.b2_mc_add_device(mc) == 0
        oks = _all_gather_obj(comm, ok)      # every device must be added before binding
        if all(oks):
            ok = lib.b2_mc_bind(mc, self.seg) == 0
            oks = _all_gather_obj(comm, ok)
        if not all(oks):
            if mc:
                lib.b2_mc_destroy(mc)
            if comm.rank == 0:
                sys.stderr.write(f"mpi4jax_b200: NVLS multicast unavailable ({native.last_error()}); "
                                 "using P2P paths only\n")
            return
        self.mc = mc
        dist.barrier(group=comm._group)

    def destroy(self) -> None:
        lib = _lib()
        if self.mc:
            lib.b2_mc_destroy(self.mc)
            self.mc = None
        if self.seg:
            lib.b2_seg_destroy(self.seg)
            self.seg = None


class NativeComm:
    """GPU side of a communicator (created collectively on first CUDA op)."""

    def __init__(self, comm: Comm):
        lib = _lib()
        setup_cuda_mpi()
        if comm.device.type != "cuda":
            raise MPIError("this process has no CUDA device; cannot communicate CUDA tensors")
        self.comm = comm
        self.device = comm.device.index
        torch.cuda.set_device(self.device)
        if lib.b2_init(self.device) != 0:
            raise MPIError(f"native init failed: {native.last_error()}")
        mode = os.environ.get("MPI4JAX_B200_HEAP", "vmm").lower()
        if mode == "vmm" and not lib.b2_vmm_supported(self.device):
            mode = "ipc"
        modes = _all_gather_obj(comm, mode)
        self.mode = "ipc" if "ipc" in modes else "vmm"
        self.want_mc = (
            self.mode == "vmm"
            and env_flag("MPI4JAX_B200_NVLS", True)
            and bool(lib.b2_multicast_supported(self.device))
            and comm.size > 1
        )
        self.want_mc = all(_all_gather_obj(comm, self.want_mc))
        devs = _all_gather_obj(comm, (socket.gethostname(), self.device))
        if len({h for h, _ in devs}) != 1:
            raise MPIError("the GPU transport needs all ranks of a communicator on one NVLink node")
        self.shared_gpu = len(set(devs)) != len(devs)   # several ranks on one GPU (testing only)
        # p2p ring slot: 16 MiB stripes give 625 GB/s on a 256 MiB sendrecv, 4 MiB ones 380 GB/s (one
        # header + credit round per 64 KiB lane stripe: profiles/r2_sweep_n8.log vs r2_p2p_n2.log).  The ring
        # area is P x 8 slots per rank -- 1 GiB at 8 ranks, 0.6 % of a B200's HBM
        slot = env_int("MPI4JAX_B200_P2P_SLOT_BYTES", 16 << 20)
        ll_cap = env_int("MPI4JAX_B200_LL_BYTES", 128 << 10)
        halo_cap = env_int("MPI4JAX_B200_HALO_BYTES", 256 << 10)
        timeout = env_float("MPI4JAX_B200_TIMEOUT", 60.0)
        ctl_bytes = int(lib.b2_layout_bytes(comm.size, slot, ll_cap, halo_cap))
        self.ctl = _Segment(comm, self.device, ctl_bytes, self.mode, want_mc=False)
        self.handle = lib.b2_comm_create(self.device, comm.rank, comm.size, self.ctl.seg,
                                         slot, ll_cap, halo_cap, timeout)
        if not self.handle:
            raise MPIError(f"native communicator creation failed: {native.last_error()}")
        # transport thresholds for THIS world size on THIS GPU model (measured table, optionally overridden by
        # a tuning file: _src/tuning.py); every rank must end up with the same numbers -- the transport
        # choice is made independently on each rank from sizes and thresholds only
        from .. import tuning

        try:
            gpu_name = torch.cuda.get_device_name(self.device)
        except Exception:                       # pragma: no cover - a name is only needed to find a table
            gpu_name = None
        self.tuning = tuning.thresholds(comm.size, gpu_name)
        seen = _all_gather_obj(comm, sorted(self.tuning.items()))
        if any(t != seen[0] for t in seen):
            raise MPIError(f"the ranks disagree on the transport thresholds (MPI4JAX_B200_TUNING_FILE?): {seen}")
        if any(self.tuning[k] != tuning.NATIVE_DEFAULTS[k] for k in ("ll_max", "oneshot_max", "nvls_min")):
            lib.b2_comm_set_tuning(self.handle, self.tuning["ll_max"], self.tuning["oneshot_max"],
                                   self.tuning["nvls_min"], 0)
        if self.tuning["bcast_mc_min"] != tuning.NATIVE_DEFAULTS["bcast_mc_min"]:
            lib.b2_comm_set_option(self.handle, b"bcast_mc_min", self.tuning["bcast_mc_min"])
        self.stage: Optional[_Segment] = None
        self._stage_half = 0
        self._retired: list = []
        self._status_pool: list = []
        self._symmetric: list = []        # (base pointer, bytes, _Segment) of symmetric_empty allocations
        self._grow_stage(_MIN_STAGE)
        if comm.size > 1:
            dist.barrier(group=comm._group)

    # -- staging ---------------------------------------------------------------
    def _grow_stage(self, total_bytes: int) -> None:
        lib = _lib()
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError(
                "mpi4jax_b200: a collective needs a larger staging buffer than is allocated, "
                "which is impossible during CUDA-graph capture. Run the function once eagerly "
                "first (mpi4jax_b200.jit does) or call mpi4jax_b200.comm_reserve(nbytes, comm=comm)."
            )
        size = _MIN_STAGE
        while size < total_bytes:
            size *= 2
        torch.cuda.synchronize()
        new = _Segment(self.comm, self.device, size, self.mode, want_mc=self.want_mc)
        lib.b2_comm_set_stage(self.handle, new.seg, new.mc)
        self._stage_half = int(lib.b2_comm_stage_half(self.handle))
        if _POISON:
            # debug mode: staging never written by a peer reads back as NaN / 0xFF.. instead of
            # stale-but-plausible data (SURVEY 5.2); the barrier keeps peers from writing early
            ptr = int(lib.b2_seg_ptr(new.seg, self.comm.rank))
            torch.as_tensor(_RawDeviceBytes(ptr, new.bytes), device=f"cuda:{self.device}").fill_(0xFF)
            torch.cuda.synchronize()
            if self.comm.size > 1:
                dist.barrier(group=self.comm._group)
        old, self.stage = self.stage, new
        if old is not None:
            # Kernels get the staging pointers BY VALUE, so a CUDA graph captured earlier keeps the old
            # segment's addresses baked into its nodes (mpi4jax_b200.jit replays them for as long as the
            # function object lives).  Unmapping here would leave them dangling on every rank; the old
            # segment therefore stays mapped until the communicator is destroyed -- the growth is
            # geometric, so the retired segments together are smaller than the live one.
            self._retired.append(old)

    def ensure_stage(self, opcode: int, blk_bytes: int) -> None:
        # same formula as b2_stage_need() (csrc/b2_collectives.cu), evaluated without leaving Python
        stride = (blk_bytes + 15) & ~15
        mult = self.comm.size if opcode in (codes.OPC_ALLTOALL, codes.OPC_SCATTER, codes.OPC_REDUCE_SCATTER) else 1
        need = stride * mult + 4096
        if need > self._stage_half:
            self._grow_stage(2 * need + 8192)

    def reserve(self, nbytes: int) -> None:
        """Make sure collectives of up to ``nbytes`` per rank (alltoall / scatter / reduce_scatter: per
        peer block times size) never have to grow the staging segment again.  Collective."""
        stride = (int(nbytes) + 15) & ~15
        need = stride * self.comm.size + 4096
        if need > self._stage_half:
            self._grow_stage(2 * need + 8192)

    @property
    def has_nvls(self) -> bool:
        return self.stage is not None and self.stage.mc is not None

    # -- plumbing ----------------------------------------------------------------
    @staticmethod
    def _stream() -> int:
        return torch.cuda.current_stream().cuda_stream

    def _check(self, rc: int, opname: str) -> None:
        if rc == 0:
            return
        msg = native.last_error()
        abort_or_raise(
            f"r{self.comm.rank} | MPI_{opname} returned error code {rc}: {msg} - aborting", rc)

    def check_device_error(self) -> None:
        buf = ctypes.create_string_buffer(512)
        code = _lib().b2_comm_check_error(self.handle, buf, 512)
        if code != 0:
            abort_or_raise(buf.value.decode(), code)

    def flush(self) -> None:
        try:
            torch.cuda.synchronize(self.device)
        except RuntimeError as exc:
            self.check_device_error()
            raise MPIError(f"CUDA failure while flushing communication: {exc}") from exc
        self.check_device_error()

    def set_tuning(self, ll_max=-1, oneshot_max=-1, nvls_min=-1, max_blocks=0) -> None:
        _lib().b2_comm_set_tuning(self.handle, ll_max, oneshot_max, nvls_min, max_blocks)

    def set_option(self, key: str, value: int) -> None:
        """Runtime switches of the native communicator: ``bcast_mc_min`` (bytes), ``nvls_pipeline`` (0/1)."""
        self._check(_lib().b2_comm_set_option(self.handle, key.encode(), int(value)), "Comm_set_option")

    def get_option(self, key: str) -> int:
        """Current value of a launch parameter: ``max_blocks``, ``sm_count``, ``bcast_mc_min``, ``nvls_pipeline``."""
        value = int(_lib().b2_comm_get_option(self.handle, key.encode()))
        if value < 0:
            raise ValueError(f"unknown communicator option {key!r}")
        return value

    @property
    def max_blocks(self) -> int:
        return self.get_option("max_blocks")

    def destroy(self) -> None:
        lib = _lib()
        try:
            torch.cuda.synchronize(self.device)
        except RuntimeError:
            pass
        if self.handle:
            lib.b2_comm_destroy(self.handle)
            self.handle = None
        if self.stage is not None:
            self.stage.destroy()
            self.stage = None
        for seg in self._retired:
            seg.destroy()
        self._retired = []
        for _, _, seg in self._symmetric:
            seg.destroy()
        self._symmetric = []
        for rec in self._status_pool:
            lib.b2_status_free(rec)
        del self._status_pool[:]
        if self.ctl is not None:
            self.ctl.destroy()
            self.ctl = None

    # -- collectives -------------------------------------------------------------
    def barrier(self) -> None:
        self._check(_lib().b2_barrier(self.handle, self._stream()), "Barrier")

    def allreduce(self, x: torch.Tensor, op_code: int, algo: int = codes.ALGO_AUTO) -> torch.Tensor:
        x, dt, op_code = _prep_reduce(x, op_code)
        out = torch.empty_like(x)
        self.ensure_stage(codes.OPC_ALLREDUCE, x.numel() * x.element_size())
        rc = _lib().b2_allreduce(self.handle, x.data_ptr(), out.data_ptr(), x.numel(), dt, op_code,
                                 algo, self._stream())
        self._check(rc, "Allreduce")
        return out

    def reduce_scatter(self, x: torch.Tensor, op_code: int, algo: int = codes.ALGO_AUTO) -> torch.Tensor:
        """MPI_Reduce_scatter_block: ``x`` is ``(size, *S)``; returns op over all ranks of block ``rank``."""
        x, dt, op_code = _prep_reduce(x, op_code)
        out = torch.empty(x.shape[1:], dtype=x.dtype, device=x.device)
        blk = out.numel()
        self.ensure_stage(codes.OPC_REDUCE_SCATTER, blk * x.element_size())
        rc = _lib().b2_reduce_scatter(self.handle, x.data_ptr(), out.data_ptr(), blk, dt, op_code, algo,
                                      self._stream())
        self._check(rc, "Reduce_scatter_block")
        return out

    # -- symmetric tensors: user memory inside the symmetric heap ---------------------------------
    def symmetric_empty(self, shape, dtype: torch.dtype) -> torch.Tensor:
        """A tensor whose storage is a symmetric segment of this communicator (same size on every rank,
        mapped into every peer and bound to an NVSwitch multicast object).  Collective.  The segment
        lives as long as the communicator."""
        shape = tuple(int(d) for d in (shape if isinstance(shape, (tuple, list, torch.Size)) else (shape,)))
        itemsize = torch.empty((), dtype=dtype).element_size()
        nbytes = max(16, itemsize * int(torch.Size(shape).numel()))
        sizes = _all_gather_obj(self.comm, nbytes)
        if len(set(sizes)) != 1:
            raise MPIError(f"symmetric_empty: every rank must ask for the same size (got {sizes} bytes)")
        torch.cuda.synchronize(self.device)
        seg = _Segment(self.comm, self.device, nbytes, self.mode, want_mc=self.want_mc)
        base = int(_lib().b2_seg_ptr(seg.seg, self.comm.rank))
        self._symmetric.append((base, seg.bytes, seg))
        raw = torch.as_tensor(_RawDeviceBytes(base, seg.bytes), device=f"cuda:{self.device}")
        return raw[: itemsize * int(torch.Size(shape).numel())].view(dtype).reshape(shape)

    def _symmetric_of(self, x: torch.Tensor):
        ptr = x.data_ptr()
        for base, nbytes, seg in self._symmetric:
            if base <= ptr and ptr + x.numel() * x.element_size() <= base + nbytes:
                return seg, ptr - base
        return None, 0

    def allreduce_inplace(self, x: torch.Tensor) -> torch.Tensor:
        """SUM-allreduce of a symmetric tensor IN PLACE, reduced inside the NVSwitch: no staging copy in,
        none out (csrc/b2_collectives.cu: b2_k_allreduce_sym)."""
        if self.comm.size == 1:
            return x
        seg, off = self._symmetric_of(x)
        if seg is None or not x.is_contiguous():
            raise ValueError("allreduce_: needs a contiguous tensor (or view) from mpi4jax_b200.symmetric_empty")
        if seg.mc is None:
            raise MPIError("allreduce_: NVLS multicast is unavailable on this communicator")
        if x.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            raise TypeError("allreduce_: the in-switch reduction supports float32, bfloat16 and float16")
        if (x.numel() * x.element_size()) % 16 or off % 16:
            raise ValueError("allreduce_: the tensor must start on a 16-byte boundary and be a multiple of 16 "
                             f"bytes long (got {x.numel() * x.element_size()} bytes at offset {off})")
        dt = codes.DTYPE_CODE[x.dtype]
        mc = int(_lib().b2_mc_ptr(seg.mc)) + off
        rc = _lib().b2_allreduce_sym(self.handle, mc, x.numel(), dt, self._stream())
        self._check(rc, "Allreduce")
        return x

    def reduce(self, x: torch.Tensor, op_code: int, root: int) -> Optional[torch.Tensor]:
        x, dt, op_code = _prep_reduce(x, op_code)
        is_root = self.comm.rank == root
        out = torch.empty_like(x) if is_root else None
        self.ensure_stage(codes.OPC_REDUCE, x.numel() * x.element_size())
        rc = _lib().b2_reduce(self.handle, x.data_ptr(), out.data_ptr() if is_root else None,
                              x.numel(), dt, op_code, root, self._stream())
        self._check(rc, "Reduce")
        return out

    def scan(self, x: torch.Tensor, op_code: int) -> torch.Tensor:
        x, dt, op_code = _prep_reduce(x, op_code)
        out = torch.empty_like(x)
        self.ensure_stage(codes.OPC_SCAN, x.numel() * x.element_size())
        rc = _lib().b2_scan(self.handle, x.data_ptr(), out.data_ptr(), x.numel(), dt, op_code,
                            self._stream())
        self._check(rc, "Scan")
        return out

    def allgather(self, x: torch.Tensor) -> torch.Tensor:
        x, lay = _layout(x)
        out = torch.empty((self.comm.size, *x.shape), dtype=x.dtype, device=x.device)
        nb = x.numel() * x.element_size()
        self.ensure_stage(codes.OPC_ALLGATHER, nb)
        self._check(_lib().b2_allgather(self.handle, x.data_ptr(), out.data_ptr(), nb, _ref(lay), self._stream()),
                    "Allgather")
        return out

    def alltoall(self, x: torch.Tensor) -> torch.Tensor:
        x, lay = _layout(x, lead=True)
        out = torch.empty(x.shape, dtype=x.dtype, device=x.device)
        nb = (x.numel() // self.comm.size) * x.element_size()
        self.ensure_stage(codes.OPC_ALLTOALL, nb)
        self._check(_lib().b2_alltoall(self.handle, x.data_ptr(), out.data_ptr(), nb, _ref(lay), self._stream()),
                    "Alltoall")
        return out

    def bcast(self, x: torch.Tensor, root: int) -> torch.Tensor:
        x = _prep(x)
        nb = x.numel() * x.element_size()
        is_root = self.comm.rank == root
        out = x if is_root else torch.empty_like(x)
        self.ensure_stage(codes.OPC_BCAST, nb)
        rc = _lib().b2_bcast(self.handle, x.data_ptr() if is_root else None,
                             None if is_root else out.data_ptr(), nb, root, None, self._stream())
        self._check(rc, "Bcast")
        return out

    def gather(self, x: torch.Tensor, root: int) -> Optional[torch.Tensor]:
        x, lay = _layout(x)
        nb = x.numel() * x.element_size()
        is_root = self.comm.rank == root
        out = (torch.empty((self.comm.size, *x.shape), dtype=x.dtype, device=x.device)
               if is_root else None)
        self.ensure_stage(codes.OPC_GATHER, nb)
        rc = _lib().b2_gather(self.handle, x.data_ptr(), out.data_ptr() if is_root else None, nb,
                              root, _ref(lay), self._stream())
        self._check(rc, "Gather")
        return out

    def scatter(self, x: torch.Tensor, root: int, out_shape, dtype) -> torch.Tensor:
        is_root = self.comm.rank == root
        out = torch.empty(out_shape, dtype=dtype, device=self.comm.device)
        nb = out.numel() * out.element_size()
        src, lay = _layout(x, lead=True) if is_root else (None, None)
        self.ensure_stage(codes.OPC_SCATTER, nb)
        rc = _lib().b2_scatter(self.handle, src.data_ptr() if is_root else None, out.data_ptr(), nb,
                               root, _ref(lay), self._stream())
        self._check(rc, "Scatter")
        return out

    # -- point to point ------------------------------------------------------------
    def _status_record(self, status: Optional[Status], itemsize: int):
        if status is None:
            return None
        rec = getattr(status, "_record", None)      # one host-mapped record per Status object
        if rec is None:
            # records of collected Status objects are reused (a Status per loop iteration must not
            # leak pinned host memory); they are freed with the communicator
            rec = self._status_pool.pop() if self._status_pool else _lib().b2_status_alloc()
            if not rec:
                raise MPIError(f"allocating a status record failed: {native.last_error()}")
            status._record = rec
            pool = self._status_pool
            weakref.finalize(status, pool.append, rec)
        return rec

    def _bind_status(self, status: Optional[Status], rec, itemsize: int) -> None:
        if status is None:
            return
        if torch.cuda.is_current_stream_capturing():
            # inside a graph the record is rewritten on every replay; read it after replay
            status._bind_native(rec, _NullEvent(self.device), itemsize)
            return
        ev = torch.cuda.Event()
        ev.record()
        status._bind_native(rec, ev, itemsize)

    def send(self, x: torch.Tensor, dest: int, tag: int) -> None:
        x = _prep(x)
        rc = _lib().b2_send(self.handle, x.data_ptr(), x.numel() * x.element_size(), dest, tag,
                            self._stream())
        self._check(rc, "Send")

    def recv(self, template: torch.Tensor, source: int, tag: int,
             status: Optional[Status]) -> torch.Tensor:
        out = torch.empty(template.shape, dtype=template.dtype, device=self.comm.device)
        rec = self._status_record(status, out.element_size())
        rc = _lib().b2_recv(self.handle, out.data_ptr(), out.numel() * out.element_size(), source, tag,
                            rec, self._stream())
        self._check(rc, "Recv")
        self._bind_status(status, rec, out.element_size())
        return out

    def sendrecv(self, sendbuf: torch.Tensor, recv_template: torch.Tensor, source: int, dest: int,
                 sendtag: int, recvtag: int, status: Optional[Status]) -> torch.Tensor:
        sendbuf = _prep(sendbuf)
        out = torch.empty(recv_template.shape, dtype=recv_template.dtype, device=self.comm.device)
        rec = self._status_record(status, out.element_size())
        rc = _lib().b2_sendrecv(self.handle, sendbuf.data_ptr(),
                                sendbuf.numel() * sendbuf.element_size(), dest, sendtag,
                                out.data_ptr(), out.numel() * out.element_size(), source, recvtag,
                                rec, self._stream())
        self._check(rc, "Sendrecv")
        self._bind_status(status, rec, out.element_size())
        return out

    # -- tensor-parallel linear: tcgen05 GEMM + in-switch allreduce (csrc/b2_gemm.cu) ----------
    def gemm_allreduce(self, x: torch.Tensor, weight: torch.Tensor) -> torch.Tensor:
        """``allreduce_SUM(x @ weight.T)`` for bf16 ``x (M, K)``, ``weight (N, K)`` in ONE kernel."""
        M, K = x.shape
        N = weight.shape[0]
        out = torch.empty((M, N), dtype=torch.bfloat16, device=x.device)
        if self.comm.size > 1:
            if not self.has_nvls:
                raise MPIError("gemm_allreduce needs NVLS multicast support")
            self.ensure_stage(codes.OPC_ALLREDUCE, M * N * 2)
        rc = _lib().b2_gemm_allreduce(self.handle, x.data_ptr(), weight.data_ptr(), out.data_ptr(), M, N, K,
                                      self._stream())
        self._check(rc, "Allreduce")
        return out

    # -- fused halo exchange ---------------------------------------------------------
    def halo_exchange(self, fields, kinds, west, east, south, north, periodic_x=True,
                      at_east_wall=False, at_north_wall=False, sw=-1, se=-1, nw=-1, ne=-1) -> None:
        """Fused single-phase 8-neighbour halo exchange (csrc/b2_halo.cu).  ``fields`` are
        float32 ``(ny, nx)`` tensors with unit inner stride and a common row pitch."""
        d = native.B2HaloDesc()
        d.nfields = len(fields)
        ny, nx = fields[0].shape
        pitch = fields[0].stride(0)
        for k, (f, kind) in enumerate(zip(fields, kinds)):
            if (f.dtype != torch.float32 or tuple(f.shape) != (ny, nx) or f.stride(1) != 1
                    or f.stride(0) != pitch):
                raise ValueError("halo_exchange needs float32 fields of one shape and row pitch")
            d.field[k] = f.data_ptr()
            d.kind[k] = {"h": 0, "u": 1, "v": 2}[kind]
        d.ny, d.nx, d.pitch = ny, nx, pitch
        d.west, d.east, d.south, d.north = west, east, south, north
        d.sw, d.se, d.nw, d.ne = sw, se, nw, ne
        d.periodic_x = int(periodic_x)
        d.at_east_wall = int(at_east_wall)
        d.at_north_wall = int(at_north_wall)
        self._check(_lib().b2_halo_exchange(self.handle, ctypes.byref(d), self._stream()), "Halo")


def _nvtx_wrap(name: str, fn):
    @functools.wraps(fn)
    def wrapped(self, *args, **kwargs):
        torch.cuda.nvtx.range_push(f"mpi4jax_b200.{name}")
        try:
            return fn(self, *args, **kwargs)
        finally:
            torch.cuda.nvtx.range_pop()

    return wrapped


#: ``MPI4JAX_B200_NVTX=1``: one NVTX range per op (visible in Nsight Systems timelines); the
#: methods are left untouched otherwise, so the fast path pays nothing (SURVEY 5.1)
NVTX_OPS = ("barrier", "allreduce", "reduce", "scan", "allgather", "alltoall", "bcast", "gather", "scatter",
            "reduce_scatter", "send", "recv", "sendrecv", "gemm_allreduce", "halo_exchange")
if env_flag("MPI4JAX_B200_NVTX", False):
    for _name in NVTX_OPS:
        setattr(NativeComm, _name, _nvtx_wrap(_name, getattr(NativeComm, _name)))


class _NullEvent:
    def __init__(self, device):
        self.device = device

    def synchronize(self):
        torch.cuda.synchronize(self.device)


def _layout(x: torch.Tensor, lead: bool = False):
    """(tensor to pass, B2Strided or None).  A non-contiguous input of a data-movement collective is
    NOT materialised by a separate torch copy kernel: its strides travel to the native kernel, which
    gathers the elements while it stages them (the fused pack of SURVEY C5).  ``lead``: dimension 0
    indexes the per-peer blocks (alltoall, scatter on the root).  Layouts the kernel cannot describe
    (more than 4 non-mergeable dimensions, overlapping / negative strides) fall back to a copy."""
    if x.numel() == 0 or (x.is_contiguous() and x.data_ptr() % 16 == 0):
        return x, None
    if x.is_contiguous():
        return x.clone(), None
    shape, stride = list(x.shape), list(x.stride())
    blk_stride = 0
    if lead:
        blk_stride = stride[0]
        shape, stride = shape[1:], stride[1:]
    dims = [(n, st) for n, st in zip(shape, stride) if n != 1]
    merged = []
    for n, st in dims:                       # merge dimensions that are contiguous with respect to each other
        if merged and merged[-1][1] == st * n:
            merged[-1] = (merged[-1][0] * n, st)
        else:
            merged.append((n, st))
    if not merged:
        merged = [(1, 1)]
    if len(merged) > 4 or any(st < 0 for _, st in merged) or blk_stride < 0:
        return x.contiguous(), None
    lay = native.B2Strided()
    lay.nd, lay.esize = len(merged), x.element_size()
    for d, (n, st) in enumerate(merged):
        lay.shape[d], lay.stride[d] = n, st
    lay.blk_stride = blk_stride
    return x, lay


def _ref(lay):
    return ctypes.byref(lay) if lay is not None else None


def _prep(x: torch.Tensor) -> torch.Tensor:
    if not x.is_contiguous():
        x = x.contiguous()
    if x.data_ptr() % 16 != 0 and x.numel() > 0:
        x = x.clone()
    return x


_BOOL_OP = {
    codes.SUM: codes.LOR, codes.MAX: codes.LOR, codes.LOR: codes.LOR, codes.BOR: codes.LOR,
    codes.PROD: codes.LAND, codes.MIN: codes.LAND, codes.LAND: codes.LAND, codes.BAND: codes.LAND,
    codes.LXOR: codes.LXOR, codes.BXOR: codes.LXOR,
}


def _prep_reduce(x: torch.Tensor, op_code: int):
    x = _prep(x)
    if x.dtype not in codes.DTYPE_CODE:
        raise TypeError(f"dtype {x.dtype} is not supported by mpi4jax_b200 reductions")
    dt = codes.DTYPE_CODE[x.dtype]
    if x.dtype == torch.bool:
        op_code = _BOOL_OP[op_code]
    elif x.dtype.is_complex and op_code not in (codes.SUM, codes.PROD):
        raise NotImplementedError("only SUM and PROD are defined for complex dtypes")
    elif x.dtype.is_floating_point and op_code not in (codes.SUM, codes.PROD, codes.MIN, codes.MAX):
        raise NotImplementedError("logical/bitwise reductions need an integer or bool dtype")
    return x, dt, op_code
